"""Static spatial adjacency stacks for the three skeleton layouts.

Mirrors the public surface of the reference generator
(`/root/reference/model/layers/graph.py:4-348`): ``Graph(layout)`` with
``get_all_adjacency() -> float64 [2, V, V]`` = (``connect``: identity + bones,
``part``: semantic left/right/limb pairs, zero diagonal), plus
``get_adjacency()`` / ``get_adjacency_type(type)``.

The reference builds the matrices from raw-skeleton joint ids and a
``use_joint`` re-indexing table; here the edges are stored directly in the
compact index space the model sees (0..V-1), which is the only form the hot
path ever consumes.  ``tests/test_layers.py`` checks every matrix against the
golden copies dumped from the reference (``tests/golden/adjacency.npz``).

Other skeletons (up to ``MAX_JOINTS`` joints) are added to the same table with
``register_layout``; every consumer of a layout name (``Graph``, the models'
``layout=`` argument, ``data.mirror``, ``DevicePrefetcher(mirror_layout=)``)
then accepts the new name.
"""
import numpy as np

# (i, j) with i < j, already in model joint order.
_EDGES = {
    "h36m": dict(
        joints=22,
        bones="0-1 0-8 1-2 2-3 4-5 4-8 5-6 6-7 8-9 8-10 9-10 9-12 9-17 10-11 12-13 13-14 14-15 "
              "14-16 17-18 18-19 19-20 19-21",
        parts="0-4 0-13 0-18 1-5 1-14 1-19 2-6 3-7 4-13 4-18 5-14 5-19 12-17 13-18 14-19 15-20 16-21",
    ),
    "cmu": dict(
        joints=25,
        bones="0-1 0-8 1-2 2-3 4-5 4-8 5-6 6-7 8-9 9-10 9-13 9-19 10-11 11-12 13-14 14-15 15-16 "
              "15-18 16-17 19-20 20-21 21-22 21-24 22-23",
        parts="0-2 0-3 0-4 0-5 0-14 0-15 0-20 0-21 1-3 1-4 1-5 1-7 1-15 1-20 2-6 4-6 4-7 4-15 4-20 "
              "4-21 5-7 5-14 5-21 13-15 13-16 13-17 13-18 13-19 13-20 14-19 14-20 14-21 15-20 15-21 "
              "16-18 16-22 17-18 17-23 18-24 19-21 19-22 19-23 19-24 22-24 23-24",
    ),
    "3dpw": dict(
        joints=23,
        bones="0-2 0-3 1-2 1-4 2-5 3-6 4-7 5-8 6-9 7-10 8-11 8-12 8-13 11-12 11-13 11-14 12-15 "
              "13-16 15-17 16-18 17-19 18-20 19-21 20-22",
        parts="0-1 0-13 0-15 1-13 1-15 3-4 3-17 3-18 4-17 4-18 6-7 6-19 6-20 7-19 7-20 9-10 12-13 "
              "15-16 17-18 19-20 21-22",
    ),
}


# the BatchNorm kernels hold the per-joint constants of a channel in one table of this many rows
MAX_JOINTS = 128


def _parse(spec):
    return [tuple(int(t) for t in e.split("-")) for e in spec.split()]


def _int(x, what):
    if isinstance(x, (bool, np.bool_)) or not isinstance(x, (int, np.integer)):
        raise TypeError(f"{what} must be an int, got {x!r}")
    return int(x)


def _edge_list(pairs, joints, what):
    out, seen = [], set()
    for e in pairs:
        if len(e) != 2:
            raise ValueError(f"{what}: {e!r} is not a pair of joint indices")
        i, j = _int(e[0], what), _int(e[1], what)
        if i == j:
            raise ValueError(f"{what}: self loop {i}-{j} (the identity is added by the graph itself)")
        if not 0 <= i < j < joints:
            raise ValueError(f"{what}: edge {i}-{j} must satisfy 0 <= i < j < joints = {joints}")
        if (i, j) in seen:
            raise ValueError(f"{what}: duplicate edge {i}-{j}")
        seen.add((i, j))
        out.append(f"{i}-{j}")
    return " ".join(out)


def register_layout(name, joints, bones, parts, mirror=None):
    """Add a skeleton layout under ``name``: ``joints`` joints (1 .. ``MAX_JOINTS``), the ``bones`` of the ``connect``
    adjacency and the semantic ``parts`` pairs, each a sequence of ``(i, j)`` with ``0 <= i < j < joints`` and no
    duplicates.  ``mirror`` is an optional ``(right, left)`` pair of equal-length, disjoint joint-index lists of the
    raw windows that ``data.mirror`` swaps; without it, mirroring the layout raises.  A name can be registered once
    and the built-in layouts cannot be replaced."""
    if not isinstance(name, str) or not name:
        raise ValueError(f"layout name must be a non-empty string, got {name!r}")
    if name in _EDGES:
        raise ValueError(f"layout {name!r} is already registered")
    joints = _int(joints, "joints")
    if not 1 <= joints <= MAX_JOINTS:
        raise ValueError(f"joints = {joints} outside 1 .. {MAX_JOINTS}")
    spec = dict(joints=joints, bones=_edge_list(bones, joints, "bones"), parts=_edge_list(parts, joints, "parts"))
    if mirror is not None:
        if len(mirror) != 2:
            raise ValueError("mirror must be a (right, left) pair of joint-index lists")
        right, left = ([_int(k, "mirror") for k in side] for side in mirror)
        if len(right) != len(left):
            raise ValueError(f"mirror: right has {len(right)} joints, left {len(left)}")
        if min(right + left, default=0) < 0:
            raise ValueError("mirror: negative joint index")
        if len(set(right)) != len(right) or len(set(left)) != len(left) or set(right) & set(left):
            raise ValueError("mirror: right and left must be disjoint lists of distinct joints")
        spec["mirror"] = (right, left)
    _EDGES[name] = spec


def mirror_lists(layout):
    """``(right, left)`` lists given to ``register_layout`` for ``layout``, or None if it was registered without."""
    return _EDGES[layout].get("mirror")


class Graph:
    """Skeleton graph of one dataset layout (``h36m`` 22 joints, ``cmu`` 25, ``3dpw`` 23, or a registered one)."""

    def __init__(self, layout="h36m"):
        if layout not in _EDGES:
            # same error class as the reference (graph.py:296-297)
            raise NotImplementedError()
        spec = _EDGES[layout]
        self.layout = layout
        self.num_joint = spec["joints"]
        self.bone_pair = [list(e) for e in _parse(spec["bones"])]
        self.part_pair = [list(e) for e in _parse(spec["parts"])]

    def _sym(self, pairs, diag):
        adj = np.eye(self.num_joint) if diag else np.zeros((self.num_joint, self.num_joint))
        for i, j in pairs:
            adj[i, j] = adj[j, i] = 1
        return adj

    def get_adjacency(self):
        return self._sym(self.bone_pair + self.part_pair, True)

    def get_adjacency_type(self, type="self"):
        if type == "self":
            return np.eye(self.num_joint)
        if type == "connect":
            return self._sym(self.bone_pair, True)
        if type == "part":
            return self._sym(self.part_pair, False)
        if type == "all":
            return self.get_adjacency()
        raise ValueError(f"Invalid graph type {type}")

    def get_all_adjacency(self):
        return np.stack([self.get_adjacency_type("connect"), self.get_adjacency_type("part")], axis=0)
