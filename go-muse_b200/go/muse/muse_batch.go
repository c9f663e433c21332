package muse

/*
#include "muse_b200.h"
*/
import "C"

import (
	"fmt"
	"runtime"
	"unsafe"
)

// Batch runs a z-normalized cross correlation between a reference series and every series of a
// comparison Group on the GPU while tracking the resulting scores (go-muse muse_batch.go:13-130).
type Batch struct {
	n           int
	ref         []float64
	batch       *C.muse_batch
	gen         uint64 // generation of the Group's device store the C batch was created on
	err         error  // what the last Run could not do (Run itself returns nil, as go-muse's does)
	Comparison  *Group
	Results     *Results
	Concurrency int
}

// Err returns the error of the last Run, or nil.  go-muse's Run cannot fail and always returns nil
// (muse_batch.go:99-130); this one can -- a CUDA error, a grouping the device store cannot key (more than 64 key
// bits) -- and keeps the signature, so a failed Run is told apart from an empty result here.
func (b *Batch) Err() error { return b.err }

// NewBatch creates a new instance with a reference timeseries, a comparison group and results.
// Errors: a comparison series of another length (muse_batch.go:24-28); a constant reference,
// "Invalid input query, Standard deviation of zero" (muse_batch.go:38-41).
func NewBatch(ref *Series, comp *Group, results *Results, cc int) (*Batch, error) {
	for _, s := range comp.series {
		if ref.Length() != s.Length() {
			return nil, fmt.Errorf("%s from comparison group series does not have the same length as the reference", s.UID())
		}
	}
	if cc < 1 {
		cc = 1
	}
	b := &Batch{ref: append([]float64(nil), ref.Values()...), Comparison: comp, Results: results, Concurrency: cc}
	// installed before anything can create the C batch: a Batch on a group that is empty now binds lazily in Run
	runtime.SetFinalizer(b, func(b *Batch) {
		if b.batch != nil {
			C.muse_batch_destroy(b.batch)
		}
	})
	if len(comp.series) == 0 {
		return b, nil
	}
	if err := b.bind(); err != nil {
		return nil, err
	}
	return b, nil
}

func (b *Batch) bind() error {
	if err := b.Comparison.syncDevice(); err != nil {
		return err
	}
	if b.batch != nil && b.gen == b.Comparison.gen {
		return nil
	}
	if b.batch != nil {
		C.muse_batch_destroy(b.batch)
		b.batch = nil
	}
	c, err := deviceContext()
	if err != nil {
		return err
	}
	rc := C.muse_batch_create(c, b.Comparison.store, (*C.double)(unsafe.Pointer(&b.ref[0])), C.int64_t(len(b.ref)), &b.batch)
	if rc != C.MUSE_OK {
		if rc == C.MUSE_ERR_STDDEV_ZERO {
			return fmt.Errorf("Invalid input query, %v", "Standard deviation of zero")
		}
		return lastError(rc)
	}
	b.gen = b.Comparison.gen
	b.n = int(C.muse_batch_fft_len(b.batch))
	return nil
}

// Run calculates the top N graphs with the highest scores; one score per distinct combination of
// the groupByLabels values, or per series when none are given.  Always returns nil, like go-muse; Err() tells
// whether the run could be carried out.
func (b *Batch) Run(groupByLabels []string) error {
	b.err = nil
	if len(b.Comparison.series) == 0 {
		return nil
	}
	if err := b.bind(); err != nil {
		b.err = err
		return nil
	}
	b.err = b.run(groupByLabels, nil, nil)
	return nil
}

// RunWhere is Run over the series of Comparison.FilterByLabelValues(labels) only, on the resident device store (no second
// store, no upload): Results end up as NewBatch(ref, <a Group of those series>, ...).Run(groupByLabels) leaves them.  When
// nothing can match -- empty labels, a key or a value no series of the group has -- it returns at once and Results are
// untouched.  Always returns nil, like Run; Err() tells whether the run could be carried out.
func (b *Batch) RunWhere(labels *Labels, groupByLabels []string) error {
	b.err = nil
	if len(b.Comparison.series) == 0 || labels == nil || labels.Len() == 0 {
		return nil
	}
	if err := b.bind(); err != nil { // uploads series added since the last call: the dictionary then knows every value
		b.err = err
		return nil
	}
	cols, ids, ok := b.Comparison.whereCols(labels)
	if !ok {
		return nil
	}
	b.err = b.run(groupByLabels, cols, ids)
	return nil
}

// run scores the bound store (whereCols / whereIDs: only the series with those label ids, muse_batch_run_where) and pushes
// the device's records through Results.Update.
func (b *Batch) run(groupByLabels []string, whereCols, whereIDs []int32) error {
	comp := b.Comparison
	r := b.Results
	cols := comp.keyCols(groupByLabels)
	topN := r.TopN
	if topN < 1 {
		return nil
	}
	scores := make([]float64, topN)
	lags := make([]int64, topN)
	idx := make([]int64, topN)
	var nOut C.int64_t
	var colPtr *C.int32_t
	if len(cols) > 0 {
		colPtr = (*C.int32_t)(unsafe.Pointer(&cols[0]))
	}
	var rc C.int
	if len(whereCols) > 0 {
		rc = C.muse_batch_run_where(b.batch, (*C.int32_t)(unsafe.Pointer(&whereCols[0])), (*C.int32_t)(unsafe.Pointer(&whereIDs[0])),
			C.int32_t(len(whereCols)), colPtr, C.int32_t(len(cols)), C.int64_t(r.MaxLag), C.int64_t(topN),
			C.double(r.Threshold), C.int32_t(r.SignFilter), C.MUSE_MODE_AUTO, 0,
			(*C.double)(unsafe.Pointer(&scores[0])), (*C.int64_t)(unsafe.Pointer(&lags[0])),
			(*C.int64_t)(unsafe.Pointer(&idx[0])), &nOut)
	} else {
		rc = C.muse_batch_run(b.batch, colPtr, C.int32_t(len(cols)), C.int64_t(r.MaxLag), C.int64_t(topN),
			C.double(r.Threshold), C.int32_t(r.SignFilter),
			(*C.double)(unsafe.Pointer(&scores[0])), (*C.int64_t)(unsafe.Pointer(&lags[0])),
			(*C.int64_t)(unsafe.Pointer(&idx[0])), &nOut)
	}
	if rc != C.MUSE_OK {
		return lastError(rc)
	}
	// the device applied the Results filter and kept the TopN best; pushing those through
	// Results.Update leaves the heap exactly as pushing every group score would
	for i := 0; i < int(nOut); i++ {
		r.Update(Score{Labels: comp.series[idx[i]].Labels(), Lag: int(lags[i]), PercentScore: scores[i]})
	}
	return nil
}
