"""Scripted episodes (ddls_b200/workload.py) in the layout the CPU oracle's batch driver takes: per episode and env-step a
template id and its mount scalars."""
import numpy as np

MOUNT_FIELDS = ('max_acceptable_jct', 'part_op_mem', 'part_dep_size', 'flow_size', 'n_mounted_workers', 'n_mounted_channels')


def script_of(wl):
    """Workload -> (template ids [B, L] int32, mount scalars [B, L] oracle MOUNT_DTYPE)."""
    from oracle.oracle import MOUNT_DTYPE
    tid = np.ascontiguousarray(wl.actions['template_id'].T, dtype=np.int32)
    mount = np.zeros(tid.shape, dtype=MOUNT_DTYPE)
    for f in MOUNT_FIELDS:
        mount[f] = wl.actions[f].T
    return tid, mount


def engine_actions(engine, tid, mount, tmap=None):
    """[B, L] script -> one ACTION_DTYPE row array per env-step; ``tmap`` maps script ids to engine template ids."""
    B, L = tid.shape
    out = []
    for s in range(L):
        a = np.zeros(B, dtype=engine.ACTION_DTYPE)
        t = tid[:, s]
        a['template_id'] = t if tmap is None else np.where(t >= 0, np.asarray(tmap, dtype=np.int32)[np.maximum(t, 0)], -1)
        for f in MOUNT_FIELDS:
            a[f] = mount[f][:, s]
        out.append(a)
    return out
