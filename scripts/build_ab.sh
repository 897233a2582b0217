#!/bin/bash
# Builds HEAD's library as madrona_b200/libmadrona_b200_A.so (git-ignored) next to
# the working tree's libmadrona_b200.so, for scripts/ab_bench.sh.
set -e
cd "$(dirname "$0")/.."
git stash -q
make -C madrona_b200 -j8 > /dev/null
cp madrona_b200/libmadrona_b200.so madrona_b200/libmadrona_b200_A.so
git stash pop -q
make -C madrona_b200 -j8 > /dev/null
ls -la madrona_b200/*.so
