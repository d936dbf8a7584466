"""Per-phase timeline of the persistent chain kernel (TT_CHAIN_TRACE=1): for every task phase, when its first task
started and its last task ended (us from the kernel's first task), the mean / max task duration, and where a task's
time goes: the mean gap before each traced event (epilogue thread 0's view; events in the order they occur).  Runs the
chain alone (pooled rows already in the workspace) and inside a whole step (pooled gather -> chain), `reps` traced
launches of each; times are means over all tasks of all launches, phase bounds medians over the launches.
GPU box only:  python scripts/chain_timeline.py [B] [P] [precision] [table] [reps]"""
import os
import subprocess
import sys

import numpy as np
import torch

os.environ["TT_CHAIN_TRACE"] = "1"
os.environ["TT_CHAIN"] = "1"
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from two_towers_overlords_b200 import TwoTowersModel, _native as N  # noqa: E402
from two_towers_overlords_b200.training import FusedTrainer  # noqa: E402

B = int(sys.argv[1]) if len(sys.argv) > 1 else 2048
P = int(sys.argv[2]) if len(sys.argv) > 2 else 512
prec = sys.argv[3] if len(sys.argv) > 3 else "bf16x3"
table = len(sys.argv) > 4 and sys.argv[4] == "table"
reps = int(sys.argv[5]) if len(sys.argv) > 5 else 5
H, Lq, Ld = 384, 32, 256
N_CTAS, SLOTS = 160, 128  # kTraceCtas, kTraceSlots (tt_step_ws.cuh)
# event kinds of tt_chain_sm100.cu (EV_*)
EVENTS = ["start", "end", "acc", "stats_in", "y_out", "y_in", "part_out", "stats_loaded", "stored", "all_in"]
NAMES = ["S", "T", "F1", "F2L", "DZ", "DX", "DW2", "DW1", "G"]

torch.manual_seed(0)
m = TwoTowersModel(projection_dim=P, precision=prec, train_table=table).cuda()
tr = FusedTrainer(m, 0.3, 1e-3, B, Lq, Ld, precision=prec, use_graph=False, ids_dtype=torch.int32,
                  mask_dtype=torch.uint8)
g = torch.Generator().manual_seed(1)
for t in tr.tok:
    if t.dtype == torch.uint8:
        t.fill_(1)
    else:
        t.copy_(torch.randint(999, 30522, t.shape, generator=g).to(t.dtype))
so = tr.step_obj
RTB, NC, NCH, NCF = (B + 127) // 128, (P + 127) // 128, (H + 127) // 128, P // 64
sms = torch.cuda.get_device_properties(0).multi_processor_count
kbt = [(B + 63) // 64, (2 * B + 63) // 64]
kcb = 8
while sum((k + kcb - 1) // kcb for k in kbt) > 48:
    kcb += 8
nch = sum((k + kcb - 1) // kcb for k in kbt)
counts = [sms, 0, 3 * RTB * NC, 3 * RTB * NCF, 3 * RTB * NC, 3 * RTB * NCH if table else 0, nch * NC * NC,
          nch * NC * NCH, sms]
offs = np.concatenate([[0], np.cumsum(counts)])


def traced(phases):
    """One traced launch -> {task: {event: us from the kernel's first event}}."""
    so.internal("trace", N_CTAS * SLOTS, 2, dtype=torch.int64).zero_()
    tr._fwd_bwd(0, phases, 0)
    torch.cuda.synchronize()
    raw = so.internal("trace", N_CTAS * SLOTS, 2, dtype=torch.int64).cpu().numpy().reshape(N_CTAS, SLOTS, 2)
    t0 = raw[:, :, 1][raw[:, :, 1] > 0].min()
    ev = {}
    for c in range(N_CTAS):
        for s in range(SLOTS):
            tag, t = int(raw[c, s, 0]), int(raw[c, s, 1])
            if t == 0:
                continue
            ev.setdefault(tag >> 4, {})[EVENTS[tag & 15]] = (t - t0) / 1e3
    return ev


def gaps(rows):
    """Mean gap before each event (from the previous event of the same task), events ordered by mean time."""
    kinds = [k for k in EVENTS if k != "start" and all(k in r for r in rows)]
    kinds.sort(key=lambda k: np.mean([r[k] - r["start"] for r in rows]))
    out, prev = [], ["start"] * len(rows)
    for k in kinds:
        d = [r[k] - r[p] for r, p in zip(rows, prev)]
        out.append(f"{k} +{np.mean(d):.1f}")
        prev = [k] * len(rows)
    return " | ".join(out)


def report(title, phases):
    for _ in range(3):
        tr._fwd_bwd(0, phases, 0)
    torch.cuda.synchronize()
    runs = [traced(phases) for _ in range(reps)]
    span = [max(r["end"] for r in ev.values() if "end" in r) for ev in runs]
    print(f"{title}: B={B} P={P} {prec} table={table}: {offs[-1]} tasks on {sms} CTAs, kcb={kcb}; {reps} traced launches, "
          f"first task start -> last task end {np.median(span):.1f} us (median; min {min(span):.1f}, max {max(span):.1f})")
    for k, nm in enumerate(NAMES):
        per_run = [[ev[i] for i in range(offs[k], offs[k + 1]) if i in ev and "start" in ev[i] and "end" in ev[i]]
                   for ev in runs]
        rows = [r for rr in per_run for r in rr]
        if not rows:
            continue
        med = lambda f: np.median([f(rr) for rr in per_run])  # noqa: E731
        dur = np.array([r["end"] - r["start"] for r in rows])
        print(f"  {nm:4s} {len(rows) // reps:4d} tasks: first start {med(lambda rr: min(r['start'] for r in rr)):6.1f}  "
              f"last start {med(lambda rr: max(r['start'] for r in rr)):6.1f}  "
              f"first end {med(lambda rr: min(r['end'] for r in rr)):6.1f}  "
              f"last end {med(lambda rr: max(r['end'] for r in rr)):6.1f}  task us mean {dur.mean():5.1f} max {dur.max():5.1f}")
        if nm == "F2L":  # the q task of a (row tile, column tile) and its p / n siblings do different work
            for role, segs in (("q", (0,)), ("p|n", (1, 2))):
                sub = [ev[i] for ev in runs for i in range(offs[k], offs[k + 1])
                       if (i - offs[k]) % 3 in segs and i in ev and "start" in ev[i] and "end" in ev[i]]
                print(f"       {role:4s} {gaps(sub)}")
        elif len(rows[0]) > 2:
            print(f"       {gaps(rows)}")


try:
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                         capture_output=True, text=True, timeout=30).stdout.strip()
except Exception:  # noqa: BLE001
    smi = torch.cuda.get_device_name(0)
print(f"device: {smi}")
tr._fwd_bwd(0, 1, 0)  # the pooled rows of slot 0, for the chain-alone launches
torch.cuda.synchronize()
report("chain alone", 2)
report("whole step (pooled gather -> chain)", 0)
