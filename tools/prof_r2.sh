# final ncu captures of the tensor-core kernels (one chunk of windows per launch), written to the directory given as $1
out=${1:?usage: tools/prof_r2.sh OUT_DIR}
mkdir -p "$out"
set -x
ncu --set full --clock-control none --import-source on -k regex:"conv_tc_kernel|cqt_ts_kernel|lognorm_split" --launch-skip 5 -c 5 -o "$out/r2_final_tc" -f python tools/profile_forward.py --reps 2 > "$out/pf.log" 2>&1
ls -la "$out" | tail -5
