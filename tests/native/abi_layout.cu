// Prints size and offset of every field of the records the kernels share with their host, and the constants they are
// built with, one line each. Built against include/simlod_abi.h by default; built with -DREFERENCE_HEADERS against the
// original project's HostDeviceInterface.h / structures.cuh it printed tests/golden/reference_abi_layout.txt, which
// tests/test_abi_and_library.py compares our output with line by line. Plain host code: nothing runs on a device.
#include <cstddef>
#include <cstdint>
#include <cstdio>
#ifdef REFERENCE_HEADERS
#include "HostDeviceInterface.h"
#include "helper_math.h"
#include "structures.cuh"
typedef Point Point_; typedef Chunk Chunk_; typedef OccupancyGrid OccupancyGrid_; typedef Node Node_;
typedef Uniforms Uniforms_; typedef Stats Stats_; typedef mat4 mat4_;
static const unsigned long long CONSTANTS[] = {MAX_POINTS_PER_NODE, POINTS_PER_CHUNK, MAX_DEPTH, GRID_NUM_CELLS / 32u, BATCH_STREAM_SIZE};
#else
#include "simlod_abi.h"
typedef SimlodPoint Point_; typedef SimlodChunk Chunk_; typedef SimlodOccupancyGrid OccupancyGrid_; typedef SimlodNode Node_;
typedef SimlodUniforms Uniforms_; typedef SimlodStats Stats_; typedef SimlodMat4 mat4_;
static const unsigned long long CONSTANTS[] = {SIMLOD_MAX_POINTS_PER_NODE, SIMLOD_POINTS_PER_CHUNK, SIMLOD_MAX_DEPTH, SIMLOD_GRID_WORDS,
                                               SIMLOD_BATCH_STREAM_SIZE};
#endif

#define SIZE(T) printf("sizeof %s %zu\n", #T, sizeof(T))
#define FIELD(T, f) printf("%s.%s %zu %zu\n", #T, #f, offsetof(T, f), sizeof(((T*)nullptr)->f))

int main() {
    const char* names[] = {"MAX_POINTS_PER_NODE", "POINTS_PER_CHUNK", "MAX_DEPTH", "GRID_WORDS", "BATCH_STREAM_SIZE"};
    for (int i = 0; i < 5; i++) printf("constant %s %llu\n", names[i], CONSTANTS[i]);
    SIZE(Point_); SIZE(Chunk_); SIZE(OccupancyGrid_); SIZE(Node_); SIZE(Uniforms_); SIZE(Stats_); SIZE(mat4_);
    FIELD(Point_, x); FIELD(Point_, y); FIELD(Point_, z); FIELD(Point_, color);
    FIELD(Chunk_, points); FIELD(Chunk_, size); FIELD(Chunk_, next);
    FIELD(OccupancyGrid_, values);
    FIELD(Node_, children); FIELD(Node_, counter); FIELD(Node_, numPoints); FIELD(Node_, level); FIELD(Node_, X); FIELD(Node_, Y);
    FIELD(Node_, Z); FIELD(Node_, countIteration); FIELD(Node_, countFlag); FIELD(Node_, name); FIELD(Node_, visible);
    FIELD(Node_, isFiltered); FIELD(Node_, isLeaf); FIELD(Node_, isLarge); FIELD(Node_, grid); FIELD(Node_, points);
    FIELD(Node_, voxelChunks); FIELD(Node_, numVoxels); FIELD(Node_, numVoxelsStored);
    FIELD(Uniforms_, width); FIELD(Uniforms_, height); FIELD(Uniforms_, time); FIELD(Uniforms_, fovy_rad); FIELD(Uniforms_, world);
    FIELD(Uniforms_, view); FIELD(Uniforms_, proj); FIELD(Uniforms_, transform); FIELD(Uniforms_, transform_updateBound);
    FIELD(Uniforms_, transformInv_updateBound); FIELD(Uniforms_, persistentBufferCapacity); FIELD(Uniforms_, momentaryBufferCapacity);
    FIELD(Uniforms_, frameCounter); FIELD(Uniforms_, boxMin); FIELD(Uniforms_, boxMax); FIELD(Uniforms_, showBoundingBox);
    FIELD(Uniforms_, showPoints); FIELD(Uniforms_, colorByNode); FIELD(Uniforms_, colorByLOD); FIELD(Uniforms_, colorWhite);
    FIELD(Uniforms_, doUpdateVisibility); FIELD(Uniforms_, doProgressive); FIELD(Uniforms_, LOD); FIELD(Uniforms_, useHighQualityShading);
    FIELD(Uniforms_, minNodeSize); FIELD(Uniforms_, pointSize); FIELD(Uniforms_, updateStats); FIELD(Uniforms_, enableEDL);
    FIELD(Uniforms_, edlStrength);
    FIELD(Stats_, frameID); FIELD(Stats_, numNodes); FIELD(Stats_, numInner); FIELD(Stats_, numLeaves); FIELD(Stats_, numNonemptyLeaves);
    FIELD(Stats_, numPoints); FIELD(Stats_, numVoxels); FIELD(Stats_, allocatedBytes_momentary); FIELD(Stats_, allocatedBytes_persistent);
    FIELD(Stats_, numVisibleNodes); FIELD(Stats_, numVisibleInner); FIELD(Stats_, numVisibleLeaves); FIELD(Stats_, numVisiblePoints);
    FIELD(Stats_, numVisibleVoxels); FIELD(Stats_, numChunksPoints); FIELD(Stats_, numChunksVoxels); FIELD(Stats_, batchletIndex);
    FIELD(Stats_, numPointsProcessed); FIELD(Stats_, numAllocatedChunks); FIELD(Stats_, chunkPoolSize); FIELD(Stats_, dbg);
    FIELD(Stats_, memCapacityReached);
    return 0;
}
