package muse

// Host-side value types of the facade: label sets, series handles, scores and the top-N collector.
// Nothing in this file touches the device.  The exported names and their behaviour are go-muse's
// (labels.go, series.go, scores.go, results.go of github.com/aouyang1/go-muse) because callers
// compile against them; the implementation is this repository's own: label sets are kept as a
// sorted pair list, the collector is a small sorted slice instead of a container/heap.

import (
	"math"
	"sort"
	"strings"
	"sync"

	"github.com/google/uuid"
)

// DefaultLabel names the label a Series receives when it is created without any.
const DefaultLabel = "uid"

// LabelMap maps label keys to label values.
type LabelMap map[string]string

type labelPair struct{ key, val string }

// Labels is an immutable label set.  Pairs are held sorted by key, so Keys() and ID() never sort
// the set itself.
type Labels struct {
	pairs []labelPair
	names []string
}

// NewLabels snapshots the map (later changes to it do not reach the set).
func NewLabels(m LabelMap) *Labels {
	ls := &Labels{pairs: make([]labelPair, 0, len(m)), names: make([]string, 0, len(m))}
	for k, v := range m {
		ls.pairs = append(ls.pairs, labelPair{k, v})
	}
	sort.Slice(ls.pairs, func(a, b int) bool { return ls.pairs[a].key < ls.pairs[b].key })
	for _, p := range ls.pairs {
		ls.names = append(ls.names, p.key)
	}
	return ls
}

// Len is the number of labels in the set.
func (ls *Labels) Len() int { return len(ls.pairs) }

// Keys lists the label keys in ascending order.  The slice is shared: do not modify it.
func (ls *Labels) Keys() []string { return ls.names }

// Get looks one key up by binary search.
func (ls *Labels) Get(key string) (string, bool) {
	i := sort.Search(len(ls.pairs), func(i int) bool { return ls.pairs[i].key >= key })
	if i < len(ls.pairs) && ls.pairs[i].key == key {
		return ls.pairs[i].val, true
	}
	return "", false
}

// ID renders "k1:v1,k2:v2" for the requested keys in ascending key order; keys the set does not
// have are skipped, no keys at all means every key.  As in go-muse the CALLER'S slice is sorted in
// place (Group.indexLabelValues relies on seeing it sorted afterwards).
func (ls Labels) ID(keys []string) string {
	if len(keys) == 0 {
		keys = ls.names
	} else if !sort.StringsAreSorted(keys) {
		sort.Strings(keys)
	}
	var sb strings.Builder
	for _, k := range keys {
		v, ok := ls.Get(k)
		if !ok {
			continue
		}
		if sb.Len() > 0 {
			sb.WriteByte(',')
		}
		sb.WriteString(k)
		sb.WriteByte(':')
		sb.WriteString(v)
	}
	return sb.String()
}

// Series is one timeseries and its label set.  The values are referenced, not copied, until the
// owning Group uploads them to the device.
type Series struct {
	vals []float64
	lab  *Labels
	uid  string
}

// NewSeries wraps y.  A nil or empty label set is replaced by {DefaultLabel: <random uuid>}.
func NewSeries(y []float64, labels *Labels) *Series {
	if labels == nil || labels.Len() == 0 {
		labels = NewLabels(LabelMap{DefaultLabel: uuid.New().String()})
	}
	return &Series{vals: y, lab: labels, uid: labels.ID(nil)}
}

// Length is the number of samples.
func (s *Series) Length() int { return len(s.vals) }

// Values exposes the samples; the facade never writes to them (Group.Roll replaces them by a new slice).
func (s *Series) Values() []float64 { return s.vals }

// Labels returns the label set given at construction.
func (s *Series) Labels() *Labels { return s.lab }

// UID identifies the series inside a Group: the ID over all of its labels.
func (s *Series) UID() string { return s.uid }

// Score is one result row; the JSON names are go-muse's wire format.
type Score struct {
	Labels       *Labels `json:"labels"`
	Lag          int     `json:"lag"`
	PercentScore float64 `json:"percentScore"`
}

func (s Score) magnitude() float64 { return math.Abs(s.PercentScore) }

// Scores is a list of Score.  The five methods below keep it usable with container/heap as a
// min-heap on |PercentScore|, which is how go-muse's callers may already hold it.
type Scores []Score

func (sc Scores) Len() int           { return len(sc) }
func (sc Scores) Less(a, b int) bool { return sc[a].magnitude() < sc[b].magnitude() }
func (sc Scores) Swap(a, b int)      { sc[a], sc[b] = sc[b], sc[a] }
func (sc *Scores) Push(v interface{}) {
	*sc = append(*sc, v.(Score))
}
func (sc *Scores) Pop() interface{} {
	last := len(*sc) - 1
	v := (*sc)[last]
	*sc = (*sc)[:last]
	return v
}

// SignFilter restricts results by the sign of the score.
type SignFilter int

// Untyped, as in go-muse, so that existing callers may also hold them in plain ints.
const (
	SignFilter_ANY = 0
	SignFilter_POS = 1
	SignFilter_NEG = -1
)

// Results collects the TopN scores by |PercentScore| among those with |Lag| <= MaxLag,
// |PercentScore| >= Threshold and the requested sign.  Safe for concurrent Update calls.  It is
// not reset between runs; Fetch empties it.
type Results struct {
	MaxLag     int
	TopN       int
	Threshold  float64
	SignFilter SignFilter

	mu   sync.Mutex
	kept Scores // ascending by magnitude; among equals the later arrival sits first
}

// NewResults builds an empty collector.
func NewResults(maxLag int, topN int, threshold float64, signFilter SignFilter) *Results {
	capHint := topN
	if capHint < 0 {
		capHint = 0
	}
	return &Results{MaxLag: maxLag, TopN: topN, Threshold: threshold, SignFilter: signFilter, kept: make(Scores, 0, capHint)}
}

func (r *Results) admits(s Score) bool {
	lag := s.Lag
	if lag < 0 {
		lag = -lag
	}
	if lag > r.MaxLag || !(s.magnitude() >= r.Threshold) { // a NaN score admits nothing
		return false
	}
	switch r.SignFilter {
	case SignFilter_ANY:
		return true
	case SignFilter_POS:
		return s.PercentScore > 0
	case SignFilter_NEG:
		return s.PercentScore < 0
	}
	return false
}

// Update offers one score.  Scores without labels are ignored.  Once TopN scores are held, a new
// one gets in only by being STRICTLY larger in magnitude than the smallest held.
func (r *Results) Update(s Score) {
	if s.Labels == nil {
		return
	}
	r.mu.Lock()
	defer r.mu.Unlock()
	if !r.admits(s) {
		return
	}
	m := s.magnitude()
	if len(r.kept) >= r.TopN {
		if r.TopN <= 0 || !(m > r.kept[0].magnitude()) {
			return
		}
		r.kept = r.kept[1:]
	}
	// first position whose magnitude is >= m: equal magnitudes already held stay behind the newcomer
	at := sort.Search(len(r.kept), func(i int) bool { return r.kept[i].magnitude() >= m })
	r.kept = append(r.kept, Score{})
	copy(r.kept[at+1:], r.kept[at:])
	r.kept[at] = s
}

// Fetch returns what is held in DESCENDING magnitude together with the mean magnitude (NaN when
// nothing is held) and leaves the collector empty.
func (r *Results) Fetch() (Scores, float64) {
	r.mu.Lock()
	defer r.mu.Unlock()
	n := len(r.kept)
	out := make(Scores, n)
	total := 0.0
	for i, s := range r.kept {
		out[n-1-i] = s
		total += s.magnitude()
	}
	r.kept = r.kept[:0]
	return out, total / float64(n)
}
