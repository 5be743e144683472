#!/bin/bash
# Burgers (main_Burgers1d.py problem) at N_domain = 16 000, N_boundary = 600 (M = 64 600), NB = 512, 8 GN steps:
# the unsharded one-GPU class path (--single) and the sharded path on 1, 2, 4, 8 GPUs (as many as the box has).
# Per-phase times are CUDA events, max over ranks (tools/dist_solve.py); GPP_TRACE adds the split of the sharded inverse
# into U = L^-T and the Theta^-1 sub-blocks, and the per-step split of the GN steps (stderr, *.trace).
# Afterwards: final loss and sol_sampled_pts of every sharded run against the one-GPU run (and the largest relative
# difference over the whole loss history, with the iteration where it occurs).
#   usage: tools/runs/r03_burgers_N16k.sh OUTDIR
set -u
OUT=${1:?output directory}
mkdir -p "$OUT"
nvidia-smi --query-gpu=index,name,power.limit,clocks.max.sm,memory.total --format=csv > "$OUT/gpus.csv"
NG=$(nvidia-smi -L | wc -l)
ARGS="--pde burgers --N 16000 --Nb 600 --NB 512 --gn_steps 8 --reps 1"
echo "GPP_TRACE=1 python tools/dist_solve.py $ARGS --single --dump-outputs $OUT/single" > "$OUT/commands.txt"
GPP_TRACE=1 python tools/dist_solve.py $ARGS --single --dump-outputs "$OUT/single" > "$OUT/single.jsonl" 2> "$OUT/single.trace"
for P in 1 2 4 8; do
  [ "$P" -le "$NG" ] || break
  CMD="python -m torch.distributed.run --nnodes=1 --nproc-per-node=$P --master-addr 127.0.0.1 --master-port 29631 tools/dist_solve.py $ARGS --dump-outputs $OUT/p$P"
  echo "GPP_TRACE=1 $CMD" >> "$OUT/commands.txt"
  GPP_TRACE=1 $CMD > "$OUT/p$P.jsonl" 2> "$OUT/p$P.trace"
done
python - "$OUT" <<'EOF'
import glob, json, os, sys
import numpy as np
out, N = sys.argv[1], 16000
band = max(1e-8, 10 * np.finfo(float).eps / 1e-5)
ref_loss = np.load(os.path.join(out, "single", "loss_hist.npy"))
ref_sol = np.load(os.path.join(out, "single", "sol.npy"))[:N]
for d in sorted(glob.glob(os.path.join(out, "p*/"))):
    loss, sol = np.load(os.path.join(d, "loss_hist.npy")), np.load(os.path.join(d, "sol.npy"))[:N]
    rel = np.abs(loss - ref_loss) / np.abs(ref_loss)
    r = dict(run=os.path.basename(d.rstrip("/")), final_loss=float(loss[-1]), final_loss_single=float(ref_loss[-1]),
             final_loss_rel=float(rel[-1]), sol_sampled_pts_rel=float(np.max(np.abs(sol - ref_sol)) / np.max(np.abs(ref_sol))),
             band=band, loss_hist_rel_max=float(rel.max()), loss_hist_rel_max_at_iter=int(rel.argmax()))
    r["final_loss_and_sol_within_band"] = r["final_loss_rel"] <= band and r["sol_sampled_pts_rel"] <= band
    print(json.dumps(r))
EOF
