package muse

/*
#include "muse_b200.h"
*/
import "C"

import (
	"fmt"
	"unsafe"
)

// RunMany scores several reference series against one comparison Group in a single call: what a loop
// of NewBatch(ref_q, comp, results_q, cc).Run(groupByLabels) computes in go-muse (muse_batch.go:23-130),
// with the store read once for up to 256 references at a time (muse_multi_run: the bounds of all of them as one
// bf16 contraction on the tensor cores).  results[q] receives the
// scores of refs[q]; a constant reference gets NewBatch's error in errs[q] and leaves results[q] untouched.
// Not part of go-muse's API: the reference builds one Batch per query.
func RunMany(refs []*Series, comp *Group, results []*Results, groupByLabels []string) (errs []error, err error) {
	return runMany(refs, comp, results, false, nil, groupByLabels)
}

// RunManyWhere is RunMany over the series of comp.FilterByLabelValues(labels) only, on the resident device store (one
// selection for every reference, no second store): results[q] ends up as RunMany on a Group of those series leaves it --
// what a loop of NewBatch(ref_q, comp, results_q, cc).RunWhere(labels, groupByLabels) computes (muse_multi_run_where).
// It makes the checks of RunMany.  When nothing can match -- empty labels, a key or a value no series of the group has --
// there is no device call: every results[q] is untouched and every errs[q] nil, as Batch.RunWhere does.
// Not part of go-muse's API.
func RunManyWhere(refs []*Series, comp *Group, results []*Results, labels *Labels, groupByLabels []string) (errs []error, err error) {
	return runMany(refs, comp, results, true, labels, groupByLabels)
}

// runMany is RunMany, or RunManyWhere when filter is set.
func runMany(refs []*Series, comp *Group, results []*Results, filter bool, labels *Labels, groupByLabels []string) (errs []error, err error) {
	if len(refs) != len(results) {
		return nil, fmt.Errorf("%d references but %d results", len(refs), len(results))
	}
	errs = make([]error, len(refs))
	if len(refs) == 0 || len(comp.series) == 0 {
		return errs, nil
	}
	n := comp.Length()
	r0 := results[0]
	rows := make([]float64, 0, len(refs)*n)
	for q, ref := range refs {
		if ref.Length() != n {
			return nil, fmt.Errorf("%s does not have the same length as the comparison group", ref.UID())
		}
		if rq := results[q]; rq.MaxLag != r0.MaxLag || rq.TopN != r0.TopN || rq.Threshold != r0.Threshold || rq.SignFilter != r0.SignFilter {
			return nil, fmt.Errorf("RunMany needs the same MaxLag, TopN, Threshold and SignFilter on every Results")
		}
		rows = append(rows, ref.Values()...)
	}
	if r0.TopN < 1 || (filter && (labels == nil || labels.Len() == 0)) {
		return errs, nil
	}
	if err := comp.syncDevice(); err != nil { // uploads series added since the last call: the dictionary then knows every value
		return nil, err
	}
	var whereCols, whereIDs []int32
	if filter {
		var ok bool
		if whereCols, whereIDs, ok = comp.whereCols(labels); !ok {
			return errs, nil
		}
	}
	c, err := deviceContext()
	if err != nil {
		return nil, err
	}
	cols := comp.keyCols(groupByLabels)
	var colPtr *C.int32_t
	if len(cols) > 0 {
		colPtr = (*C.int32_t)(unsafe.Pointer(&cols[0]))
	}
	topN := r0.TopN
	scores := make([]float64, len(refs)*topN)
	lags := make([]int64, len(refs)*topN)
	idx := make([]int64, len(refs)*topN)
	nOut := make([]int64, len(refs))
	var rc C.int
	if filter {
		rc = C.muse_multi_run_where(c, comp.store, (*C.double)(unsafe.Pointer(&rows[0])), C.int64_t(len(refs)), C.int64_t(n),
			(*C.int32_t)(unsafe.Pointer(&whereCols[0])), (*C.int32_t)(unsafe.Pointer(&whereIDs[0])), C.int32_t(len(whereCols)),
			colPtr, C.int32_t(len(cols)), C.int64_t(r0.MaxLag), C.int64_t(topN), C.double(r0.Threshold),
			C.int32_t(r0.SignFilter), C.MUSE_MODE_AUTO,
			(*C.double)(unsafe.Pointer(&scores[0])), (*C.int64_t)(unsafe.Pointer(&lags[0])),
			(*C.int64_t)(unsafe.Pointer(&idx[0])), (*C.int64_t)(unsafe.Pointer(&nOut[0])))
	} else {
		rc = C.muse_multi_run(c, comp.store, (*C.double)(unsafe.Pointer(&rows[0])), C.int64_t(len(refs)), C.int64_t(n),
			colPtr, C.int32_t(len(cols)), C.int64_t(r0.MaxLag), C.int64_t(topN), C.double(r0.Threshold),
			C.int32_t(r0.SignFilter), C.MUSE_MODE_AUTO,
			(*C.double)(unsafe.Pointer(&scores[0])), (*C.int64_t)(unsafe.Pointer(&lags[0])),
			(*C.int64_t)(unsafe.Pointer(&idx[0])), (*C.int64_t)(unsafe.Pointer(&nOut[0])))
	}
	if rc != C.MUSE_OK {
		return nil, lastError(rc)
	}
	for q := range refs {
		if nOut[q] < 0 {
			errs[q] = fmt.Errorf("Invalid input query, %v", "Standard deviation of zero")
			continue
		}
		for i := 0; i < int(nOut[q]); i++ {
			k := q*topN + i
			results[q].Update(Score{Labels: comp.series[idx[k]].Labels(), Lag: int(lags[k]), PercentScore: scores[k]})
		}
	}
	return errs, nil
}
