#!/bin/sh
# Link-compatibility check ("existing callers link unchanged"): compile the reference's OWN tutorial
# tutorials/minimal/minimal.cpp, untouched and against the reference's OWN headers, and link it against
# libembree4_b200.so instead of libembree4.so.  Only the resulting binaries are kept, in oracle/_ref/link_compat with the
# other reference build products (git-ignored); no reference source enters the repo.  Runs only where the reference exists;
# elsewhere the binaries built before are used (tests/test_link_compat.py).  Our host drivers are in tests/link_compat/.
set -e
cd "$(dirname "$0")"
REF=${EMBREE_REFERENCE:-/root/reference}
GEN=_ref/gen_rel/include/embree4
[ -f "$REF/tutorials/minimal/minimal.cpp" ] && [ -d "$GEN" ] || { echo "reference not present: keeping prebuilt binary"; exit 0; }
# -lembree4 resolves to libembree4_b200.so through this alias; the binaries record the library's soname
# (libembree4_b200.so) and find it through their rpath, $ORIGIN/../../../embree_b200/csrc
OUT=_ref/link_compat
HOST=../tests/link_compat
GOLD=../tests/golden
mkdir -p $OUT
ln -sf ../../../embree_b200/csrc/libembree4_b200.so $OUT/libembree4.so
g++ -O1 -std=c++11 -I"$REF/include" -I"$GEN" -o $OUT/embree_minimal "$REF/tutorials/minimal/minimal.cpp" \
    -L$OUT -lembree4 -Wl,-rpath,'$ORIGIN/../../../embree_b200/csrc'
echo built oracle/_ref/link_compat/embree_minimal

# BASELINE configs[0]: the reference's tutorial device code tutorials/triangle_geometry/triangle_geometry_device.cpp (cube +
# ground plane, rtcTraversableIntersect1 + rtcTraversableOccluded1 per pixel in its own tile loop), compiled untouched
# together with the reference's sys / tasking sources it needs and OUR small host driver (tutorial_host.cpp: what
# tutorial.cpp would provide), linked (a) against libembree4_b200.so -> oracle/_ref/link_compat/embree_triangle_geometry (runs on the GPU
# box) and (b) against the unmodified reference library -> the golden frame tests/golden/triangle_geometry_160x120.raw.
GENR=_ref/gen_rel
INC="-I$REF -I$REF/include -I$GENR/include -I$GENR/include/embree4 -I$GENR -DTASKING_INTERNAL"
SYS="$REF/common/sys/sysinfo.cpp $REF/common/sys/alloc.cpp $REF/common/sys/thread.cpp $REF/common/sys/mutex.cpp $REF/common/sys/condition.cpp
     $REF/common/sys/barrier.cpp $REF/common/sys/estring.cpp $REF/common/sys/regression.cpp $REF/common/tasking/taskschedulerinternal.cpp
     $REF/common/math/constants.cpp $REF/tutorials/common/alloc/alloc.cpp"
if [ ! -x $OUT/embree_triangle_geometry ] || [ $HOST/tutorial_host.cpp -nt $OUT/embree_triangle_geometry ]; then
  g++ -O1 -std=c++17 -w $INC -o $OUT/embree_triangle_geometry $HOST/tutorial_host.cpp "$REF/tutorials/triangle_geometry/triangle_geometry_device.cpp" $SYS \
      -L$OUT -lembree4 -lpthread -Wl,-rpath,'$ORIGIN/../../../embree_b200/csrc'
  echo built oracle/_ref/link_compat/embree_triangle_geometry
fi
if [ -f _ref/libembree4.so.4 ] && [ ! -f $GOLD/triangle_geometry_160x120.raw ]; then
  g++ -O1 -std=c++17 -w $INC -o $OUT/ref_triangle_geometry $HOST/tutorial_host.cpp "$REF/tutorials/triangle_geometry/triangle_geometry_device.cpp" $SYS \
      -L_ref -l:libembree4.so.4 -lpthread -Wl,-rpath,'$ORIGIN/..'
  $OUT/ref_triangle_geometry $GOLD/triangle_geometry_160x120.raw 160 120 4
  rm -f $OUT/ref_triangle_geometry
fi

# BASELINE configs[3]a: the reference's tutorial device code tutorials/hair_geometry/hair_geometry_device.cpp (hair sets converted with
# rtcSetGeometryTessellationRate / rtcSetGeometryEnableFilterFunctionFromArguments, per pixel a path of rtcTraversableIntersect1 and
# rtcTraversableOccluded1 with its transparency-accumulating occlusion filter), compiled untouched with OUR host driver hair_host.cpp
# (procedural fur ball: round linear / flat Bezier / round Bezier hair), linked (a) against libembree4_b200.so ->
# oracle/_ref/link_compat/embree_hair_geometry and (b) against the unmodified reference -> golden frames tests/golden/hair_geometry_<type>_96x72.raw.
if [ ! -x $OUT/embree_hair_geometry ] || [ $HOST/hair_host.cpp -nt $OUT/embree_hair_geometry ]; then
  g++ -O1 -std=c++17 -w $INC -o $OUT/embree_hair_geometry $HOST/hair_host.cpp "$REF/tutorials/hair_geometry/hair_geometry_device.cpp" $SYS \
      -L$OUT -lembree4 -lpthread -Wl,-rpath,'$ORIGIN/../../../embree_b200/csrc'
  echo built oracle/_ref/link_compat/embree_hair_geometry
fi
if [ -f _ref/libembree4.so.4 ] && [ ! -f $GOLD/hair_geometry_2_96x72.raw ]; then
  g++ -O1 -std=c++17 -w $INC -o $OUT/ref_hair_geometry $HOST/hair_host.cpp "$REF/tutorials/hair_geometry/hair_geometry_device.cpp" $SYS \
      -L_ref -l:libembree4.so.4 -lpthread -Wl,-rpath,'$ORIGIN/..'
  for t in 0 1 2; do $OUT/ref_hair_geometry $GOLD/hair_geometry_${t}_96x72.raw 96 72 4 $t 3000; done
  rm -f $OUT/ref_hair_geometry
fi

# BASELINE configs[3]b: the reference's tutorial device code tutorials/dynamic_scene/dynamic_scene_device.cpp (DYNAMIC | ROBUST scene of a plane
# and 20 spheres with per-geometry build qualities, all vertices rewritten and re-committed every frame), compiled untouched with OUR host
# driver dynamic_host.cpp, linked (a) against libembree4_b200.so -> oracle/_ref/link_compat/embree_dynamic_scene and (b) against the unmodified reference ->
# golden frames tests/golden/dynamic_scene_160x120_<frame>.raw.
if [ ! -x $OUT/embree_dynamic_scene ] || [ $HOST/dynamic_host.cpp -nt $OUT/embree_dynamic_scene ]; then
  g++ -O1 -std=c++17 -w $INC -o $OUT/embree_dynamic_scene $HOST/dynamic_host.cpp "$REF/tutorials/dynamic_scene/dynamic_scene_device.cpp" $SYS \
      -L$OUT -lembree4 -lpthread -Wl,-rpath,'$ORIGIN/../../../embree_b200/csrc'
  echo built oracle/_ref/link_compat/embree_dynamic_scene
fi
if [ -f _ref/libembree4.so.4 ] && [ ! -f $GOLD/dynamic_scene_160x120_2.raw ]; then
  g++ -O1 -std=c++17 -w $INC -o $OUT/ref_dynamic_scene $HOST/dynamic_host.cpp "$REF/tutorials/dynamic_scene/dynamic_scene_device.cpp" $SYS \
      -L_ref -l:libembree4.so.4 -lpthread -Wl,-rpath,'$ORIGIN/..'
  $OUT/ref_dynamic_scene $GOLD/dynamic_scene_160x120 160 120 4 3
  rm -f $OUT/ref_dynamic_scene
fi

# Point primitives: the reference's tutorial device code tutorials/point_geometry/point_geometry_device.cpp (three sets of 512 sphere /
# disc / oriented-disc points over a ground plane, closest hit + shadow ray per pixel), compiled untouched with tutorial_host.cpp (camera of
# point_geometry.cpp:23-24), linked (a) against libembree4_b200.so -> oracle/_ref/link_compat/embree_point_geometry and (b) against the unmodified reference ->
# the golden frame tests/golden/point_geometry_160x120.raw.
PCAM="-DCAMERA_FROM=0.0f,2.0f,7.0f"
if [ ! -x $OUT/embree_point_geometry ] || [ $HOST/tutorial_host.cpp -nt $OUT/embree_point_geometry ]; then
  g++ -O1 -std=c++17 -w $INC $PCAM -o $OUT/embree_point_geometry $HOST/tutorial_host.cpp "$REF/tutorials/point_geometry/point_geometry_device.cpp" $SYS \
      -L$OUT -lembree4 -lpthread -Wl,-rpath,'$ORIGIN/../../../embree_b200/csrc'
  echo built oracle/_ref/link_compat/embree_point_geometry
fi
if [ -f _ref/libembree4.so.4 ] && [ ! -f $GOLD/point_geometry_160x120.raw ]; then
  g++ -O1 -std=c++17 -w $INC $PCAM -o $OUT/ref_point_geometry $HOST/tutorial_host.cpp "$REF/tutorials/point_geometry/point_geometry_device.cpp" $SYS \
      -L_ref -l:libembree4.so.4 -lpthread -Wl,-rpath,'$ORIGIN/..'
  $OUT/ref_point_geometry $GOLD/point_geometry_160x120.raw 160 120 4
  rm -f $OUT/ref_point_geometry
fi
