# builds the library of the CURRENT csrc/ into variants/<name>.so (experiments: several builds timed in one GPU visit, tools/gpu_variants.sh);
# sources and flags are agarcl_b200/build.py's, $EXTRA adds nvcc flags
set -eo pipefail
cd "$(dirname "$0")/.."
mkdir -p variants
python -c 'import shlex, subprocess, sys; sys.path.insert(0, "agarcl_b200"); import build
subprocess.check_call(build.nvcc_command(sys.argv[1], shlex.split(sys.argv[2]), verbose=True))' "variants/$1.so" "${EXTRA:-}" 2>&1 \
  | grep -A2 "k_stepENS\|error" | grep "stack\|Used\|error"
