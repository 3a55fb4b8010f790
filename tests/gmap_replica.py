"""A plain-Python restatement of the GPU-resident keypoint map (csrc/gmap.cu), for tests.

It follows the oracle's Map (src/mymap.cpp, src/keypoint.cpp:23-32, updateMap) and adds what the oracle does not keep:
the update that wrote each entry (its tag), the export order and the storable-position rule.  Every float operation is a
numpy float32 operation, so it rounds as the fp32 device code does (no FMA).

- position: R p + T as ((r0 x + r1 y) + r2 z) + t, then createKeypoint's int(trunc(v / 10)) * 10;
- block: getBlockID, int(roundf(v / 10000)) * 10000 per axis (half away from zero), 21 bits each;
- admission: rejected when an entry of the block lies within 800 mm and is at least as salient (<=); otherwise an entry at
  the same lattice position is overwritten in place (it takes the new update's tag), else the keypoint is appended;
- blocks in creation order, entries of a block in insertion order;
- a position is storable when every transformed, unsnapped coordinate is finite and within +-STORABLE_MM; other
  keypoints are skipped, and they are not dropped ones.
"""
import math

import numpy as np

f32 = np.float32
PREC = 10000
LATTICE = f32(10.0)
REJECT_MM = f32(800.0)
STORABLE_MM = f32(2.1e9)


def roundf(v):
    """C roundf of a float32: half away from zero"""
    v = float(v)
    return int(math.copysign(math.floor(abs(v) + 0.5), v))


def snap(v):
    """Keypoint::createKeypoint: int(trunc(v / 10)) * 10"""
    return f32(int(math.trunc(float(f32(v) / LATTICE))) * 10)


def block_coord(v):
    return roundf(f32(v) / f32(PREC))


def block_id(x, y, z):
    key = 0
    for v in (x, y, z):
        key = (key << 21) | ((block_coord(v) * PREC) & 0x1FFFFF)
    return key


def transform(xyz, pose):
    """R p + T in fp32 with the map update's rounding; pose = row-major 3 x 4 (None = identity)"""
    xyz = np.asarray(xyz, f32).reshape(-1, 3)
    if pose is None:
        return xyz.copy()
    P = np.asarray(pose, f32).reshape(3, 4)
    x, y, z = xyz[:, 0], xyz[:, 1], xyz[:, 2]
    with np.errstate(invalid="ignore", over="ignore"):
        return np.stack([((P[r, 0] * x + P[r, 1] * y) + P[r, 2] * z) + P[r, 3] for r in range(3)], axis=1).astype(f32)


def storable(xyz):
    with np.errstate(invalid="ignore"):
        return np.all(np.abs(np.asarray(xyz, f32)) <= STORABLE_MM, axis=-1)


class Map:
    """blocks: block id -> list of entries [x, y, z, ratio, desc (6,) uint64, tag]"""

    def __init__(self):
        self.blocks = {}
        self.updates = 0

    def __len__(self):
        return sum(len(b) for b in self.blocks.values())

    def add(self, xyz, ratio, desc, pose=None):
        """one map update (bshot_gmap_add): every keypoint in order.  Returns the number of keypoints skipped as not storable"""
        w = transform(xyz, pose)
        ratio = np.asarray(ratio, f32).reshape(-1)
        desc = np.asarray(desc, np.uint64).reshape(-1, 6)
        if len(w) == 0:
            return 0
        tag, skipped = self.updates, 0
        ok = storable(w)
        for i in range(len(w)):
            if not ok[i]:
                skipped += 1
                continue
            e = [snap(w[i, 0]), snap(w[i, 1]), snap(w[i, 2]), ratio[i], desc[i].copy(), tag]
            blk = self.blocks.setdefault(block_id(e[0], e[1], e[2]), [])
            reject, same = False, None
            for k, q in enumerate(blk):
                dx, dy, dz = e[0] - q[0], e[1] - q[1], e[2] - q[2]
                if np.sqrt((dx * dx + dy * dy) + dz * dz) < REJECT_MM and e[3] <= q[3]:
                    reject = True
                if same is None and (q[0], q[1], q[2]) == (e[0], e[1], e[2]):
                    same = k
            if reject:
                continue
            if same is None:
                blk.append(e)
            else:
                blk[same] = e
        self.updates += 1
        return skipped

    def _cube(self, pos, rng):
        pos = np.asarray(pos, f32).reshape(3)
        rng = f32(rng)
        return [(roundf((pos[a] - rng) / f32(PREC)), roundf((pos[a] + rng) / f32(PREC))) for a in range(3)]

    def probes(self, pos, rng):
        """blocks getKeypoints visits around pos"""
        c = self._cube(pos, rng)
        return max(0, c[0][1] - c[0][0] + 1) * max(0, c[1][1] - c[1][0] + 1) * max(0, c[2][1] - c[2][0] + 1)

    def get(self, pos, rng):
        """Map::getKeypoints: entries of the blocks of the +-rng cube, x outermost, z innermost -> (xyz, desc, tags)"""
        (x0, x1), (y0, y1), (z0, z1) = self._cube(pos, rng)
        out = []
        for bx in range(x0, x1 + 1):
            for by in range(y0, y1 + 1):
                for bz in range(z0, z1 + 1):
                    out += self.blocks.get(block_id(f32(bx * PREC), f32(by * PREC), f32(bz * PREC)), [])
        return _arrays(out)

    def export(self):
        """gmap_export's map order: blocks in ascending lattice coordinates -> (xyzr, desc, tags)"""
        out = []
        for blk in sorted((b for b in self.blocks.values() if b), key=lambda b: tuple(block_coord(v) for v in b[0][:3])):
            out += blk
        xyz, desc, tags = _arrays(out)
        ratio = np.array([e[3] for e in out], f32).reshape(-1, 1)
        return np.concatenate([xyz, ratio], axis=1), desc, tags


def _arrays(entries):
    xyz = np.array([e[:3] for e in entries], f32).reshape(-1, 3)
    desc = np.array([e[4] for e in entries], np.uint64).reshape(-1, 6)
    tags = np.array([e[5] for e in entries], np.uint32)
    return xyz, desc, tags
