"""Reading and writing the committed fixtures of tests/golden.

A fixture stores what a computation returned, kept small:
  * inputs are not stored: they are drawn again from their seeds here (`intree_inputs`, `nll_analysis_inputs`) and
    checked against the SHA-256 the fixture recorded of the arrays the computation was given;
  * volumes the tests compare with a tolerance are stored on a fixed, seeded sample of their voxels (`Fixture.sample`
    takes the same sample of a computed volume); volumes compared bit for bit are stored whole;
  * an array identical to an earlier one is stored once.
"""
import hashlib
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
N_SAMPLE = 4096

# v1_tta.npz / v1_notta.npz: which part of the 182x218x182 result each entry holds; the argmax is stored as packed
# bits on the voxels of `v1_seg_sample`
V1_LATTICE = np.s_[::6, ::6, ::6]          # class-1 probability on a stride-6 lattice
V1_BLOCK = np.s_[68:100, 88:120, 68:100]   # both probabilities, dense 32^3 block


def digest(a) -> str:
    a = np.ascontiguousarray(a)
    return hashlib.sha256(("%s %s " % (a.dtype.str, a.shape)).encode() + a.tobytes()).hexdigest()


def v1_seg_sample(shape):
    """A seeded half of the voxels.  Planes or lattices would follow the stride-2 structure of the network's output
    (the no-TTA foreground fraction is 0.591 over the volume, 0.604 over even z planes)."""
    return np.random.default_rng(0).random(shape, dtype=np.float32) < 0.5


def save_v1(path, seg, probs, **extra):
    m = v1_seg_sample(seg.shape)
    np.savez_compressed(path, seg_bits=np.packbits(seg[m]), shape=np.array(seg.shape), seg_sample_sha256=np.array(digest(m)),
                        p1_lattice=probs[1][V1_LATTICE].astype(np.float32), p1_block=probs[1][V1_BLOCK].astype(np.float32),
                        p0_block=probs[0][V1_BLOCK].astype(np.float32), fg_frac=np.array([seg[m].mean()]), **extra)


def load_v1(path):
    """-> dict of the stored arrays plus `seg_sample` (boolean volume) and `seg` (the argmax on those voxels)."""
    g = dict(np.load(path))
    m = v1_seg_sample(tuple(int(s) for s in g["shape"]))
    assert digest(m) == str(g["seg_sample_sha256"]), "the seeded voxel sample differs from the one the fixture stores"
    g["seg_sample"], g["seg"] = m, np.unpackbits(g["seg_bits"])[: int(m.sum())]
    return g


class Fixture(dict):
    def __init__(self, arrays, index, shape):
        super().__init__(arrays)
        self._index, self._shape = index, shape

    def sample(self, a):
        """The stored voxel sample of a volume of the fixture's shape."""
        a = np.asarray(a)
        assert a.shape == self._shape, (a.shape, self._shape)
        return a.reshape(-1)[self._index]


def save(path, arrays, inputs, sampled, seed=0):
    """arrays: name -> array to store; inputs: name -> array as the computation saw it (digest only); sampled: names of
    volumes stored on the voxel sample (all of one shape)."""
    shape = {np.shape(arrays[k]) for k in sampled}
    assert len(shape) == 1, shape
    shape = shape.pop()
    index = np.sort(np.random.default_rng(seed).choice(int(np.prod(shape)), size=N_SAMPLE, replace=False)).astype(np.int32)
    out = {"sample_index": index, "sample_shape": np.array(shape),
           "input_names": np.array(sorted(inputs)), "input_sha256": np.array([digest(inputs[k]) for k in sorted(inputs)])}
    seen = {digest(v): k for k, v in inputs.items()}
    alias_names, alias_targets = [], []
    for k, v in arrays.items():
        v = np.asarray(v)
        d = digest(v)
        if v.size > 64 and d in seen and (k in sampled or seen[d] not in sampled):
            alias_names.append(k); alias_targets.append(seen[d])
            continue
        seen.setdefault(d, k)
        out[k] = v.reshape(-1)[index] if k in sampled else v
    out["alias_names"], out["alias_targets"] = np.array(alias_names, dtype=str), np.array(alias_targets, dtype=str)
    out["sampled_names"] = np.array(sorted(sampled))
    np.savez_compressed(path, **out)


def load(path, inputs) -> Fixture:
    """Stored arrays plus the regenerated inputs (each checked against its recorded digest); aliases resolved, sampled
    names already sampled."""
    f = np.load(path)
    index, shape = f["sample_index"], tuple(int(s) for s in f["sample_shape"])
    arrays = {k: f[k] for k in f.files}
    for name, d in zip(f["input_names"].tolist(), f["input_sha256"].tolist()):
        assert digest(inputs[name]) == d, "regenerated input %s differs from the one the fixture was made from" % name
        arrays[name] = inputs[name]
    sampled = set(f["sampled_names"].tolist())
    for name, target in zip(f["alias_names"].tolist(), f["alias_targets"].tolist()):
        a = arrays[target]
        arrays[name] = a.reshape(-1)[index] if name in sampled and target not in sampled else a
    return Fixture(arrays, index, shape)


def intree() -> Fixture:
    return load(os.path.join(HERE, "intree_v1.npz"), intree_inputs())


def nll_analysis() -> Fixture:
    return load(os.path.join(HERE, "nll_analysis_v1.npz"), nll_analysis_inputs())


# ------------------------------------------------------------------------------------------------
# seeded inputs
# ------------------------------------------------------------------------------------------------
def stage1_inputs(seed=7, shape=(40, 46, 38), k=5):
    """Seeded stage-1 inputs: a target, k registered references, a rough brain mask, a valid-score mask."""
    rng = np.random.default_rng(seed)
    g = np.stack(np.meshgrid(*[np.linspace(-1, 1, s) for s in shape], indexing="ij"))
    brain = ((g ** 2).sum(0) < 0.8).astype("float32")
    base = (100 + 30 * g[0] + 20 * np.sin(3 * g[1]) * g[2]).astype("float32")
    refs = [(base * rng.uniform(0.8, 1.2) + rng.normal(0, 8, shape)).astype("float32") * brain for _ in range(k)]
    target = (base + rng.normal(0, 8, shape)).astype("float32")
    target[12:16, 20:25, 15:19] += 80.0                          # a hyper-intense lesion
    target *= brain
    valid = (brain * (rng.random(shape) > 0.1)).astype("float32")
    return target, refs, brain, valid


def masked_z_score(x, mask):
    """z-score over mask > 0 with numpy.ma statistics: bit for bit what the reference's z_score returned on the
    fixture's volumes, as float32 (its digest in intree_v1.npz checks this)."""
    m = np.ma.masked_array(x, mask=1 - mask)
    return ((x - m.mean()) / max(m.std(), 0.00001)).astype(np.float32)


def intree_inputs():
    """Everything intree_v1.npz's computations were given, in the order make_golden_intree.py draws it."""
    target, refs, brain, valid = stage1_inputs()
    rng = np.random.default_rng(11)
    sparks = (rng.random((30, 34, 28)) > 0.8).astype("float32")
    shape = (33, 40, 29)
    xs = [np.clip(rng.normal(0.5, 0.35, size=shape), 0, 1).astype(np.float32) for _ in range(5)]
    xs[2][:4] = 0.5
    m = (rng.random(shape) > 0.3).astype(np.float32)
    a = (rng.random((20, 20, 20)) > 0.6).astype("float32")
    b = (rng.random((20, 20, 20)) > 0.6).astype("float32")
    rng2 = np.random.default_rng(31)
    gm = [(rng2.random(target.shape) > 0.35).astype("float32") for _ in refs]
    for x in gm:
        x[5:9] = 0                                               # a slab no reference covers -> NaN
    speck = valid.copy()
    speck[2:4, 3:6, 4:6] = 1.0                                   # sparks outside the brain, to be filtered away
    speck[36:39, 40:43, 30:34] = 1.0
    zt = masked_z_score(target, brain)
    return {"in_target": target, "in_refs": np.stack(refs), "in_brain": brain, "in_valid": valid, "sparks_in": sparks,
            "ens_x": np.stack(xs), "ens_mask": m, "dice_in": np.stack([a, b]), "gmask": np.stack(gm), "cf_in": speck,
            "z_target": zt, "zscore_masked": zt, "z_refs": np.stack([masked_z_score(r, brain) for r in refs])}


def nll_analysis_inputs():
    """The case nll_analysis_v1.npz's run was given: target, k references, their brain masks and tissue labels."""
    rng = np.random.default_rng(23)
    shape, k = (44, 52, 40), 6
    g = np.stack(np.meshgrid(*[np.linspace(-1, 1, s) for s in shape], indexing="ij"))
    r2 = (g ** 2).sum(0)
    base = (100 + 25 * g[0] + 15 * np.cos(2 * g[1]) * g[2]).astype("float32")
    brains, tissues, refs = [], [], []
    for i in range(k):
        rad = 0.78 + 0.04 * rng.random()
        brain = (r2 < rad).astype("float32")
        # tissue labels 0..3 (background / cerebrum / cerebellum + brainstem / cortex), slightly different per reference
        t = np.zeros(shape, "float32")
        t[r2 < rad] = 3
        t[r2 < rad - 0.12] = 1
        t[(r2 < rad - 0.05) & (g[2] < -0.35 + 0.03 * rng.random()) & (g[1] < 0.1)] = 2
        img = ((base * rng.uniform(0.85, 1.15) + rng.normal(0, 7, shape)) * brain).astype("float32")
        refs.append(img); brains.append(brain); tissues.append(t)
    target = (base + rng.normal(0, 7, shape)).astype("float32")
    target[14:18, 22:27, 20:24] += 70.0                              # lesion in the cerebrum
    target[20:23, 12:15, 6:9] += 60.0                                # lesion in the cerebellum (median-filtered region)
    target *= (r2 < 0.8)
    return {"in_target": target, "in_refs": np.stack(refs), "in_label1": np.stack(brains),
            "in_label2": np.stack(tissues).astype(np.uint8)}
