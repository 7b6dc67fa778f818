// bridge.go — the thin cgo layer between the reference's Go package `core` and the B200
// library (include/rs_knn.h -> librs_knn_b200.so).  This file is what a maintainer of
// Oneaccount1/recommend-sys adds; it could not be compiled in the build image (no Go
// toolchain), so every behaviour it relies on is exercised through the same C ABI by the
// Python mirror (recommend-sys_b200/core.py) and the C++ mirror (host/core.hpp).
//
// cgo rules honoured here:
//   - C never retains a Go pointer: every slice is borrowed for the duration of one call
//     (rs_knn_fit / rs_knn_predict_batch copy to the device before returning);
//   - goroutines migrate between OS threads, so the library binds the CUDA device on every
//     entry (api.cu: enter());
//   - Go `int` is 64-bit: inner ids are narrowed to int32 when marshalled;
//   - the handle lives in an UNEXPORTED field so gob (core/dump.go:11-43, used by Copy in
//     core/eval.go:29-30) neither serialises nor aliases it.
package core

/*
#cgo CFLAGS: -I${SRCDIR}/../../../include
#cgo LDFLAGS: -L${SRCDIR}/../.. -lrs_knn_b200 -Wl,-rpath,${SRCDIR}/../..
#include <stdlib.h>
#include "rs_knn.h"
*/
import "C"

import (
	"fmt"
	"reflect"
	"runtime"
	"unsafe"
)

// simEnum maps a Sim func value to the library's enum by comparing code pointers
// (core/sim.go:7 makes Sim a plain func type; the device cannot call back into Go).
// Any other function is an error: there is no CPU fallback.
func simEnum(s Sim) C.int32_t {
	p := reflect.ValueOf(s).Pointer()
	switch p {
	case reflect.ValueOf(Cosine).Pointer():
		return C.RS_SIM_COSINE
	case reflect.ValueOf(MSD).Pointer():
		return C.RS_SIM_MSD
	case reflect.ValueOf(Pearson).Pointer():
		return C.RS_SIM_PEARSON
	case reflect.ValueOf(PearsonBaseline).Pointer():
		return C.RS_SIM_PEARSON_BASELINE
	}
	panic("core: the CUDA KNN supports the built-in similarities only (Cosine, MSD, Pearson, PearsonBaseline)")
}

func knnTypeEnum(t string) C.int32_t {
	switch t {
	case basic:
		return C.RS_KNN_BASIC
	case centered:
		return C.RS_KNN_CENTERED
	case zScore:
		return C.RS_KNN_ZSCORE
	case baseline:
		return C.RS_KNN_BASELINE
	}
	panic("core: unknown KNN type " + t)
}

// check panics on a non-zero status: the reference has no error returns on this path
// (core/base.go:68-74 panics, core/base.go:26-54 type assertions panic).
func check(rc C.int32_t) {
	if rc != C.RS_OK {
		panic(fmt.Sprintf("rs_knn error %d: %s", int(rc), C.GoString(C.rs_last_error())))
	}
}

type deviceKNN struct{ h *C.rs_knn }

func newDeviceKNN(p Parameters, knnType string) *deviceKNN {
	var cp C.rs_knn_params
	check(C.rs_knn_params_default(&cp))
	cp.sim = simEnum(p.GetSim("sim", MSD))
	cp.knn_type = knnTypeEnum(knnType)
	cp.k = C.int32_t(p.GetInt("k", 40))
	cp.min_k = C.int32_t(p.GetInt("mink", 1))
	cp.device = C.int32_t(p.GetInt("device", -1))
	if p.GetString("pearsonMode", "exact") == "sums" {
		cp.pearson_mode = C.RS_PEARSON_SUMS
	}
	switch p.GetString("simPath", "auto") {
	case "tensor":
		cp.sim_path = C.RS_PATH_TENSOR
	case "stream":
		cp.sim_path = C.RS_PATH_STREAM
	}
	if p.GetString("store", "matrix") == "topk" {
		cp.store = C.RS_STORE_TOPK
	}
	cp.topk = C.int32_t(p.GetInt("topk", p.GetInt("k", 40)))
	cp.row_begin = C.int64_t(p.GetInt("rowBegin", 0))
	cp.row_end = C.int64_t(p.GetInt("rowEnd", 0))
	cp.shrinkage = C.double(p.GetFloat64("shrinkage", 0))
	// sharding over the GPUs of one box (rs_knn.h: symmetric slabs for RS_STORE_TOPK, cyclic row
	// shards for RS_STORE_MATRIX); 0 = this handle computes everything
	cp.shard_count = C.int32_t(p.GetInt("shardCount", 0))
	cp.shard_index = C.int32_t(p.GetInt("shardIndex", 0))
	d := &deviceKNN{}
	check(C.rs_knn_create(&cp, &d.h))
	runtime.SetFinalizer(d, func(d *deviceKNN) { d.close() })
	return d
}

func (d *deviceKNN) close() {
	if d.h != nil {
		C.rs_knn_destroy(d.h)
		d.h = nil
	}
}

func i32(p []int32) *C.int32_t {
	if len(p) == 0 {
		return nil
	}
	return (*C.int32_t)(unsafe.Pointer(&p[0]))
}

func f64(p []float64) *C.double {
	if len(p) == 0 {
		return nil
	}
	return (*C.double)(unsafe.Pointer(&p[0]))
}

func (d *deviceKNN) fit(left, right []int32, rating []float64, nLeft, nRight int, globalMean float64,
	leftBias, rightBias []float64, globalBias float64) {
	check(C.rs_knn_fit(d.h, i32(left), i32(right), f64(rating), C.int64_t(len(rating)),
		C.int32_t(nLeft), C.int32_t(nRight), C.double(globalMean), f64(leftBias), f64(rightBias),
		C.double(globalBias)))
	runtime.KeepAlive(left)
	runtime.KeepAlive(right)
	runtime.KeepAlive(rating)
}

// update adds ratings (inner ids, in call order) to the fitted model: it becomes the Fit of the union (rs_knn_update).
func (d *deviceKNN) update(left, right []int32, rating []float64, nLeft, nRight int, globalMean float64) {
	check(C.rs_knn_update(d.h, i32(left), i32(right), f64(rating), C.int64_t(len(rating)), C.int32_t(nLeft),
		C.int32_t(nRight), C.double(globalMean)))
	runtime.KeepAlive(left)
	runtime.KeepAlive(right)
	runtime.KeepAlive(rating)
}

// baselineALS is the EXTENSION behind Parameters["baseline"] = "als" (BASELINE.json config 3): ALS
// baseline estimates computed on the device instead of BaseLine.Fit's sequential SGD
// (core/base.go:135-163).  Returns (userBias, itemBias); the global bias is the global mean.
func baselineALS(device int, users, items []int32, rating []float64, nUsers, nItems int, globalMean,
	regU, regI float64, nEpochs int) ([]float64, []float64) {
	ub, ib := make([]float64, nUsers), make([]float64, nItems)
	check(C.rs_baseline_als(C.int32_t(device), i32(users), i32(items), f64(rating), C.int64_t(len(rating)),
		C.int32_t(nUsers), C.int32_t(nItems), C.double(globalMean), C.double(regU), C.double(regI),
		C.int32_t(nEpochs), f64(ub), f64(ib)))
	return ub, ib
}

// setK forwards Parameters["k"] / ["mink"], which the reference reads at Predict time
// (core/knn.go:80-81), to a fitted handle.
func (d *deviceKNN) setK(k, minK int) { check(C.rs_knn_set_k(d.h, C.int32_t(k), C.int32_t(minK))) }

// Cyclic row shards (one estimator per GPU, Parameters["shardCount"] >= 2 with the matrix kept):
// peerExport returns the 64-byte CUDA IPC handle + offset of this shard's matrix, peerImport
// attaches all shards' matrices (gathered by whatever transport joins the processes), mirror pulls
// the triangle this shard did not compute over NVLink.  With all shards in ONE process
// (goroutine per GPU, like the reference's nJobs) peerImportLocal takes the handles directly.
func (d *deviceKNN) peerExport() ([64]byte, int64) {
	var hb [64]byte
	var off C.int64_t
	check(C.rs_knn_peer_export(d.h, (*C.uchar)(unsafe.Pointer(&hb[0])), &off))
	return hb, int64(off)
}

func (d *deviceKNN) peerImport(handles [][64]byte, offsets []int64) {
	flat := make([]byte, 64*len(handles))
	for i := range handles {
		copy(flat[64*i:], handles[i][:])
	}
	check(C.rs_knn_peer_import(d.h, C.int32_t(len(handles)), (*C.uchar)(unsafe.Pointer(&flat[0])),
		(*C.int64_t)(unsafe.Pointer(&offsets[0]))))
}

func (d *deviceKNN) peerImportLocal(peers []*deviceKNN) {
	hs := make([]*C.rs_knn, len(peers))
	for i, p := range peers {
		hs[i] = p.h
	}
	check(C.rs_knn_peer_import_local(d.h, C.int32_t(len(hs)), &hs[0]))
}

func (d *deviceKNN) mirror() { check(C.rs_knn_mirror(d.h)) }

// predictBatchShardedDevice: every shard gets the FULL test set (device pointers), answers the pairs whose left
// row it owns and leaves +0.0 elsewhere (a cold-start pair is answered by shard index % shardCount); an int64 SUM
// all-reduce of the bit patterns over the shards (NCCL) then holds the complete prediction vector on every GPU.
func (d *deviceKNN) predictBatchShardedDevice(dLeft, dRight unsafe.Pointer, n int, dOut unsafe.Pointer) {
	check(C.rs_knn_predict_batch_sharded_device(d.h, (*C.int32_t)(dLeft), (*C.int32_t)(dRight), C.int64_t(n),
		(*C.double)(dOut)))
}

// recommendShardedDevice: every shard gets the same queries (device pointers) and writes its PARTIAL lists
// ids[n][nTop] / scores[n][nTop]: the targets it owns for right queries, the whole list of the left queries whose row
// it owns.  All-gather them and unite them with rs_knn_topk_union_device (groups of at most 2048 / nTop lists).
func (d *deviceKNN) recommendShardedDevice(side int, dQueries unsafe.Pointer, n, nTop int, dIDs, dScores unsafe.Pointer) {
	check(C.rs_knn_recommend_sharded_device(d.h, C.int32_t(side), (*C.int32_t)(dQueries), C.int64_t(n), C.int32_t(nTop),
		(*C.int32_t)(dIDs), (*C.double)(dScores)))
}

// scoreAllShardedDevice: the score rows out[n][nTargets] of this shard, +0.0 in the cells it does not answer; an
// int64 SUM all-reduce of the bit patterns over the shards assembles rs_knn_score_all.
func (d *deviceKNN) scoreAllShardedDevice(side int, dQueries unsafe.Pointer, n int, dOut unsafe.Pointer) {
	check(C.rs_knn_score_all_sharded_device(d.h, C.int32_t(side), (*C.int32_t)(dQueries), C.int64_t(n),
		(*C.double)(dOut)))
}

func (d *deviceKNN) predictBatch(left, right []int32) []float64 {
	out := make([]float64, len(left))
	check(C.rs_knn_predict_batch(d.h, i32(left), i32(right), C.int64_t(len(left)), f64(out)))
	return out
}

// Query sides of rs_knn_recommend (enum rs_side).
const (
	sideLeft  = 0
	sideRight = 1
)

// recommend: ids / scores are [len(queries)][nTop], row-major.
func (d *deviceKNN) recommend(side int, queries []int32, nTop int) ([]int32, []float64) {
	ids := make([]int32, len(queries)*nTop)
	scores := make([]float64, len(queries)*nTop)
	if len(queries) == 0 {
		return ids, scores
	}
	check(C.rs_knn_recommend(d.h, C.int32_t(side), i32(queries), C.int64_t(len(queries)), C.int32_t(nTop), i32(ids),
		f64(scores)))
	return ids, scores
}

// recommendGiven: queries given as rating lists — list b is ids[ptr[b]:ptr[b+1]] (inner ids of the target side) with
// ratings vals[...], in the caller's order (rs_knn_recommend_given).  ids / scores are [len(ptr)-1][nTop], row-major.
func (d *deviceKNN) recommendGiven(side int, ptr []int64, ids []int32, vals []float64, nTop int) ([]int32, []float64) {
	n := len(ptr) - 1
	outIDs := make([]int32, n*nTop)
	outScores := make([]float64, n*nTop)
	if n <= 0 {
		return outIDs, outScores
	}
	if len(ids) == 0 { // every list empty: the library still wants valid pointers
		ids, vals = []int32{0}, []float64{0}
	}
	check(C.rs_knn_recommend_given(d.h, C.int32_t(side), (*C.int64_t)(unsafe.Pointer(&ptr[0])), i32(ids), f64(vals),
		C.int64_t(n), C.int32_t(nTop), i32(outIDs), f64(outScores)))
	return outIDs, outScores
}

// pinnedInt32 / pinnedFloat64: page-locked host memory of the library's per-process cache (rs_knn_host_alloc) viewed
// as a Go slice, for callers that stage large batches themselves: copies from and to such memory run at full PCIe
// speed.  The memory is C memory (no Go pointers in it); release returns the block to the cache.
func pinnedInt32(n int) (s []int32, release func()) {
	var p unsafe.Pointer
	check(C.rs_knn_host_alloc(C.size_t(n*4), &p))
	return unsafe.Slice((*int32)(p), n), func() { C.rs_knn_host_free(p) }
}

func pinnedFloat64(n int) (s []float64, release func()) {
	var p unsafe.Pointer
	check(C.rs_knn_host_alloc(C.size_t(n*8), &p))
	return unsafe.Slice((*float64)(p), n), func() { C.rs_knn_host_free(p) }
}

func (d *deviceKNN) simsRows(row0, nrows, n int) []float64 {
	out := make([]float64, nrows*n)
	check(C.rs_knn_sims_rows(d.h, C.int64_t(row0), C.int64_t(nrows), f64(out)))
	return out
}

func (d *deviceKNN) topK(k, rows int) ([]int32, []float64) {
	idx := make([]int32, rows*k)
	sim := make([]float64, rows*k)
	check(C.rs_knn_topk(d.h, C.int32_t(k), i32(idx), f64(sim)))
	return idx, sim
}

func (d *deviceKNN) means(n int) []float64 {
	out := make([]float64, n)
	check(C.rs_knn_means(d.h, f64(out)))
	return out
}

func (d *deviceKNN) stddevs(n int) []float64 {
	out := make([]float64, n)
	check(C.rs_knn_stddevs(d.h, f64(out)))
	return out
}
