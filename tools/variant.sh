# Build a variant of one translation unit with extra -D flags into libmcmcn_<name>.so (same ABI; A/B with tools/ab.sh):
#   bash tools/variant.sh <name> -DMCMCN_DEBUG_BOUNDS                     (the tcgen05 step kernel, mcmcn_sets_tc.cu)
#   UNIT=mcmcn_sets_logit bash tools/variant.sh <name> -DMY_SWITCH=1 ...   (a switch added to the source for the A/B)
set -e
name=$1; shift
unit=${UNIT:-mcmcn_sets_tc}
root=$(cd "$(dirname "$0")/.." && pwd)
csrc=$root/mcmc-for-nested-data_b200/csrc
/usr/local/cuda/bin/nvcc -gencode arch=compute_100a,code=sm_100a -lineinfo -O3 -std=c++17 -I $root/include -I $csrc -Xcompiler -fPIC "$@" \
  -c $csrc/$unit.cu -o /tmp/${unit}_$name.o
objs=$(ls $csrc/build/*.o | grep -v $unit.o)
/usr/local/cuda/bin/nvcc -shared --cudart shared -o $root/mcmc-for-nested-data_b200/libmcmcn_$name.so $objs /tmp/${unit}_$name.o -ldl
echo built libmcmcn_$name.so
