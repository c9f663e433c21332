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

// Sharded comparison groups: one process per GPU of a box (MUSE_DEVICE = local rank), each holding a contiguous
// block of the group's series; the reference is given to every process.  go-muse has no such mode -- its Batch.Run
// walks one in-memory Group (muse_batch.go:99-130) -- so this file is an addition, not a mirror: the scores,
// the group max before the filter (muse_batch.go:87-89), the filter (results.go:46-52) and the top-N
// (results.go:54-87) of the WHOLE group come out of every process identical to a single-process Run.
//
// A step is one call, Batch.RunSharded: the kernels that produce a shard's records store them into every process's
// receive buffer over NVLink peer memory and the merge runs on the device (muse_batch_run_exchange_ex); there is no
// collective library underneath.  Setup needs one out-of-band exchange of 64 bytes per process (Handle /
// OpenPeers), e.g. over the launcher's rendezvous.

// ExchangeHandleBytes is the size of the handle every process publishes to its peers.
const ExchangeHandleBytes = 64

// Exchange is this process's end of the peer-memory exchange.
type Exchange struct {
	x     *C.muse_exchange
	rank  int
	world int
}

// NewExchange creates the receive buffers for `capacity` records per peer and step: at least TopN for runs without
// groupByLabels, at least the number of label groups a shard can hold for grouped runs.
func NewExchange(rank, world, capacity int) (*Exchange, error) {
	c, err := deviceContext()
	if err != nil {
		return nil, err
	}
	if world < 1 || rank < 0 || rank >= world {
		return nil, fmt.Errorf("muse_b200: rank %d of %d", rank, world)
	}
	e := &Exchange{rank: rank, world: world}
	if rc := C.muse_exchange_create(c, C.int32_t(rank), C.int32_t(world), C.int64_t(capacity), &e.x); rc != C.MUSE_OK {
		return nil, lastError(rc)
	}
	runtime.SetFinalizer(e, func(e *Exchange) { e.Close() })
	return e, nil
}

// Handle returns the 64 bytes the other processes need to map this process's receive buffers.
func (e *Exchange) Handle() ([]byte, error) {
	h := make([]byte, ExchangeHandleBytes)
	if rc := C.muse_exchange_ipc_handle(e.x, unsafe.Pointer(&h[0])); rc != C.MUSE_OK {
		return nil, lastError(rc)
	}
	return h, nil
}

// OpenPeers maps every process's buffers; handles[r] is what rank r's Handle returned.
func (e *Exchange) OpenPeers(handles [][]byte) error {
	if len(handles) != e.world {
		return fmt.Errorf("muse_b200: %d handles for %d ranks", len(handles), e.world)
	}
	all := make([]byte, 0, e.world*ExchangeHandleBytes)
	for r, h := range handles {
		if len(h) != ExchangeHandleBytes {
			return fmt.Errorf("muse_b200: handle of rank %d has %d bytes", r, len(h))
		}
		all = append(all, h...)
	}
	if rc := C.muse_exchange_open_peers(e.x, unsafe.Pointer(&all[0])); rc != C.MUSE_OK {
		return lastError(rc)
	}
	return nil
}

// Close releases the buffers (peers must have stopped stepping).
func (e *Exchange) Close() {
	if e.x != nil {
		C.muse_exchange_destroy(e.x)
		e.x = nil
	}
}

// SetShard declares this Group to be the block of a sharded group that starts at series index `first` of the whole,
// and fixes the label dictionary: for every label key the complete list of its values, IDENTICAL on every
// process, so that the int32 ids the device groups by mean the same labels everywhere.  Call before the first
// NewBatch on the group.
func (g *Group) SetShard(first int64, dictionary map[string][]string) {
	g.sharded = true
	g.shardFirst = first
	g.fixedDict = dictionary
	if g.store != nil { // re-encode with the fixed ids
		C.muse_group_destroy(g.store)
		g.store = nil
		g.uploaded = 0
	}
}

// ShardScore is one score of the whole sharded group.  Index counts series over all shards in rank order; Labels is
// set when that series lives in this process's shard (the other processes hold the rest).
type ShardScore struct {
	Index        int64
	Lag          int
	PercentScore float64
	Labels       *Labels
}

// RunSharded is Batch.Run over the whole sharded group: every process calls it the same number of times with the same
// groupByLabels and Results settings, and every process gets the same scores back, best first (results.go:54-87).
func (b *Batch) RunSharded(e *Exchange, groupByLabels []string) ([]ShardScore, error) {
	comp := b.Comparison
	if len(comp.series) == 0 {
		return nil, errNoSeries
	}
	if err := b.bind(); err != nil {
		return nil, err
	}
	r := b.Results
	if r.TopN < 1 {
		return nil, nil
	}
	cols := comp.keyCols(groupByLabels)
	scores := make([]float64, r.TopN)
	lags := make([]int64, r.TopN)
	idx := make([]int64, r.TopN)
	var nOut C.int64_t
	var colPtr *C.int32_t
	if len(cols) > 0 {
		colPtr = (*C.int32_t)(unsafe.Pointer(&cols[0]))
	}
	rc := C.muse_batch_run_exchange_ex(b.batch, e.x, colPtr, C.int32_t(len(cols)), C.int64_t(r.MaxLag), C.int64_t(r.TopN),
		C.double(r.Threshold), C.int32_t(r.SignFilter), C.MUSE_MODE_AUTO,
		(*C.double)(unsafe.Pointer(&scores[0])), (*C.int64_t)(unsafe.Pointer(&lags[0])),
		(*C.int64_t)(unsafe.Pointer(&idx[0])), &nOut)
	if rc != C.MUSE_OK {
		return nil, lastError(rc)
	}
	out := make([]ShardScore, int(nOut))
	for i := range out {
		out[i] = ShardScore{Index: idx[i], Lag: int(lags[i]), PercentScore: scores[i]}
		if local := idx[i] - comp.shardFirst; local >= 0 && local < int64(len(comp.series)) {
			out[i].Labels = comp.series[local].Labels()
		}
	}
	return out, nil
}

// RunManySharded is RunMany over the whole sharded group (without groupByLabels): refs[q] is scored against the series of
// every process, and scores[q] -- identical on every process, best first, filled as RunSharded fills its result -- is what a
// single-process RunMany over the whole group puts into results[q].  results supply the settings (the same MaxLag, TopN,
// Threshold and SignFilter on every Results) and are left untouched.  A constant reference gets NewBatch's error in errs[q].
// Every process calls it with the same references and settings; a process whose shard holds no series takes part all the
// same.  One call runs the queries in steps of up to 256, each one exchange step (muse_multi_run_exchange).
func RunManySharded(e *Exchange, refs []*Series, comp *Group, results []*Results) (errs []error, scores [][]ShardScore, err error) {
	if len(refs) != len(results) {
		return nil, nil, fmt.Errorf("%d references but %d results", len(refs), len(results))
	}
	errs = make([]error, len(refs))
	scores = make([][]ShardScore, len(refs))
	if len(refs) == 0 {
		return errs, scores, nil
	}
	if len(comp.series) == 0 && comp.n == 0 { // an empty shard: its store takes the references' length
		comp.n = refs[0].Length()
	}
	n := comp.Length()
	r0 := results[0]
	rows := make([]float64, 0, len(refs)*n)
	for q, ref := range refs {
		if ref.Length() != n {
			return nil, nil, fmt.Errorf("%s does not have the same length as the comparison group", ref.UID())
		}
		if rq := results[q]; rq.MaxLag != r0.MaxLag || rq.TopN != r0.TopN || rq.Threshold != r0.Threshold || rq.SignFilter != r0.SignFilter {
			return nil, nil, fmt.Errorf("RunManySharded needs the same MaxLag, TopN, Threshold and SignFilter on every Results")
		}
		rows = append(rows, ref.Values()...)
	}
	if r0.TopN < 1 {
		return errs, scores, nil
	}
	if err := comp.syncDevice(); err != nil {
		return nil, nil, err
	}
	topN := r0.TopN
	sc := make([]float64, len(refs)*topN)
	lags := make([]int64, len(refs)*topN)
	idx := make([]int64, len(refs)*topN)
	nOut := make([]int64, len(refs))
	rc := C.muse_multi_run_exchange(comp.store, e.x, (*C.double)(unsafe.Pointer(&rows[0])), C.int64_t(len(refs)), C.int64_t(n),
		C.int64_t(r0.MaxLag), C.int64_t(topN), C.double(r0.Threshold), C.int32_t(r0.SignFilter), C.MUSE_MODE_AUTO,
		(*C.double)(unsafe.Pointer(&sc[0])), (*C.int64_t)(unsafe.Pointer(&lags[0])),
		(*C.int64_t)(unsafe.Pointer(&idx[0])), (*C.int64_t)(unsafe.Pointer(&nOut[0])))
	if rc != C.MUSE_OK {
		return nil, nil, lastError(rc)
	}
	for q := range refs {
		if nOut[q] < 0 {
			errs[q] = fmt.Errorf("Invalid input query, %v", "Standard deviation of zero")
			continue
		}
		out := make([]ShardScore, int(nOut[q]))
		for i := range out {
			k := q*topN + i
			out[i] = ShardScore{Index: idx[k], Lag: int(lags[k]), PercentScore: sc[k]}
			if local := idx[k] - comp.shardFirst; local >= 0 && local < int64(len(comp.series)) {
				out[i].Labels = comp.series[local].Labels()
			}
		}
		scores[q] = out
	}
	return errs, scores, nil
}
